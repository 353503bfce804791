"""--no-pairing (MM_F_INDEPEND_SEG, worker_for map.c:458-498): the two reads of a pair are flipped per pe_ori as for a joint
pair, then each is mapped on its own, and the records still print as a pair.  So the exact oracle is this build's own
single-segment path: mate 1 must map as mm_map_frag(n_segs=1) of mate 1 under its own name, mate 2 as mm_map_frag(n_segs=1)
of revcomp(mate 2) with qs/qe/rev flipped back, and no hit may carry proper_frag.  The CLI's records must equal those of the
single-end runs on r1 and on revcomp(r2) once the pairing fields are set aside."""
import ctypes as C
import hashlib
import os
import subprocess
import numpy as np
import pytest
import _libs as L
from test_gpu_api import Reg1, StepHead, _hit
from test_gpu_paths import data  # noqa: F401  (fixture: repeat family, overlapping mates, z-drop cuts)

pytestmark = pytest.mark.gpu
SYN = os.path.join(L.ROOT, "build", "mmsynth")
NEW = os.path.join(L.ROOT, "build", "minimap2-b200")
MM_F_CIGAR, MM_F_OUT_SAM, MM_F_FRAG_MODE, MM_F_INDEPEND_SEG = 0x004, 0x008, 0x2000, 0x20000

# size and sha256 of the --no-pairing CLI outputs of test_cli_equals_single_end, for machines without oracle/_ref/minimap2_B
# source: this project's output on a B200, recorded where no reference build was available; the test also holds every record,
# field by field, to the single-end runs, so these guard against regressions rather than prove parity with the reference
CLI_DIGESTS = {
    "--no-pairing -ax sr -t 8 ref.fa r1.fq r2.fq":
        {"bytes": 3415672, "sha256": "e597f5bc51c8bc8ec501de0eb0390c2f0f8a91bf8f12bab4191c00e084493803"},
    "--no-pairing -ax sr --secondary=yes -t 8 ref.fa r1.fq r2.fq":
        {"bytes": 4040679, "sha256": "4c573c789dffcefb219dd066f138e3f168be933fba8f4338931dc07d1fbda962"},
    "--no-pairing -ax sr --cs --MD -t 8 ref.fa r1.fq r2.fq":
        {"bytes": 3518525, "sha256": "65c979d8ce51ef8e8dc54c2620e9c6af1536001984feb28155006f9c9bd90d7e"},
    "--no-pairing -cx sr -t 8 ref.fa r1.fq r2.fq":
        {"bytes": 1184499, "sha256": "85c5ece5959f203a869a4480b3f84c6fb22db94067480a3c6d2a5f81d221c968"},
}


def _fastq(name, seq, qual=None):
    return b"@" + name + b"\n" + seq + b"\n+\n" + (qual if qual is not None else b"I" * len(seq)) + b"\n"


def _read_fq(fn):
    ls = open(fn, "rb").read().split(b"\n")
    return [(ls[i][1:].split()[0], ls[i + 1], ls[i + 3]) for i in range(0, len(ls) - 3, 4)]


def _write_rc(src, dst):
    """the reads of src reverse-complemented (qualities reversed), names kept"""
    with open(dst, "wb") as f:
        for n, s, q in _read_fq(src):
            f.write(_fastq(n, L.revcomp(s), q[::-1]))


# ---------------------------------------------------------------------------------------------------- device layer

def test_device_flips_from_table():
    """mmg_batch_t.flip: single-read fragments whose flips come from a table chain exactly as the same reads uploaded
    already reverse-complemented (K1-K3 and the re-chain pass see one-segment units)."""
    import airlift_b200.api as api
    from test_oracle_vs_ref import _mk_ref, _frags
    rng = np.random.default_rng(11)
    refseqs = _mk_ref(rng, n_ctg=2, ln=60000)
    ctx = api.Context(0)
    idx = api.Index(ctx, refseqs, 11, 21)
    try:
        mapped = _frags(rng, refseqs, 300, True)  # [m1, revcomp(m2)]
        opt = api.sr_opt()
        units = [[s] for f in mapped for s in (f[0], L.revcomp(f[1]))]      # the reads as read, one per unit
        flips = np.array([j for _ in mapped for j in (0, 1)], dtype=np.uint8)
        want_b, keep_w = api.Context.make_batch([[s] for f in mapped for s in f])
        want = api.chains_to_py(ctx.seed_chain_batch(idx, opt, want_b))
        got_b, keep_g = api.Context.make_batch(units)
        ctx.batch_upload(opt, got_b, flips)
        got = api.chains_to_py(ctx.seed_chain_resident(idx, opt, True))
        for k in ("n_u", "n_a", "rep_len", "n_mini", "rechained", "u_off", "a_off", "mini_off"):
            assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k
        assert np.asarray(got["u"]).tobytes() == np.asarray(want["u"]).tobytes()
        assert np.asarray(got["a"]).tobytes() == np.asarray(want["a"]).tobytes()
        assert np.array_equal(got["mini_pos"], want["mini_pos"])
        assert int(np.asarray(want["n_u"]).sum()) > 300
        with pytest.raises(ValueError):
            ctx.batch_upload(opt, got_b, flips[:-1])
    finally:
        idx.close()
        ctx.close()


# ---------------------------------------------------------------------------------------------------- library API

class Api:
    def __init__(self, ref, preset):
        import bench
        self.bench = bench
        lib = self.lib = bench.load_lib()
        lib.mm_map_frag.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.c_int),
                                    C.POINTER(C.POINTER(Reg1)), C.c_void_p, C.POINTER(bench.MapOptFull), C.c_char_p]
        lib.mm_tbuf_init.restype = C.c_void_p
        lib.mm_tbuf_destroy.argtypes = [C.c_void_p]
        self.ipt, self.opt = bench.IdxOpt(), bench.MapOptFull()
        lib.mm_set_opt(None, C.byref(self.ipt), C.byref(self.opt))
        lib.mm_set_opt(preset, C.byref(self.ipt), C.byref(self.opt))
        self.opt.flag |= MM_F_CIGAR | MM_F_OUT_SAM
        rd = lib.mm_idx_reader_open(str(ref).encode(), C.byref(self.ipt), None)
        self.mi = lib.mm_idx_reader_read(rd, 4)
        lib.mm_idx_reader_close(rd)
        lib.mm_mapopt_update(C.byref(self.opt), self.mi)
        self.tb = lib.mm_tbuf_init()

    def opt_with(self, flag):
        o = self.bench.MapOptFull()
        C.memmove(C.byref(o), C.byref(self.opt), C.sizeof(o))
        o.flag |= flag
        return o

    def read_batch(self, fns, opt):
        arr = (C.c_char_p * len(fns))(*[str(f).encode() for f in fns])
        reader = self.lib.mm_b200_open_reads(len(fns), arr)
        b = self.lib.mm_b200_read_batch(reader, C.byref(opt), 10**9)
        self.lib.mm_b200_close_reads(reader)
        return b

    @staticmethod
    def batch_hits(b):
        """{read: ([hit tuple + proper_frag], rep_len)} of a mapped batch"""
        h = C.cast(b, C.POINTER(StepHead)).contents
        return [([_hit(h.reg[r][i]) + (h.reg[r][i].bits >> 13 & 1,) for i in range(h.n_reg[r])], h.rep_len[r]) for r in range(h.n_seq)]

    def map_frag(self, name, seqs, opt, flip_qlen=None):
        n = len(seqs)
        arr = (C.c_char_p * n)(*seqs)
        qlens = (C.c_int * n)(*[len(s) for s in seqs])
        n_regs = (C.c_int * n)()
        regs = (C.POINTER(Reg1) * n)()
        self.lib.mm_map_frag(self.mi, n, qlens, arr, n_regs, regs, self.tb, C.byref(opt), name)
        out = [[_hit(regs[j][i], flip_qlen) + (regs[j][i].bits >> 13 & 1,) for i in range(n_regs[j])] for j in range(n)]
        rep_len = C.cast(self.tb, C.POINTER(C.c_int))[0]  # mm_tbuf_t: {rep_len, frag_gap}
        return out, rep_len

    def close(self):
        self.lib.mm_tbuf_destroy(self.tb)
        self.lib.mm_idx_destroy(self.mi)


def _check_independent(api, r1, r2, flip2, every=1):
    """map r1/r2 as pairs with MM_F_INDEPEND_SEG through mm_b200_map_batch; every `every`-th pair must equal
    mm_map_frag(n_segs=1) of each mate (mate 2 reverse-complemented when flip2, its hits flipped back).  Returns the batch hits,
    the number of hits checked and the path counters of the batch call."""
    opt = api.opt_with(MM_F_INDEPEND_SEG)
    b = api.read_batch([r1, r2], opt)
    pc = (C.c_uint64 * 8)()
    api.lib.mm_b200_path_counts(api.mi, pc, 1)
    assert api.lib.mm_b200_map_batch(api.mi, C.byref(opt), 8, b, 0) == 0
    api.lib.mm_b200_path_counts(api.mi, pc, 1)
    got = api.batch_hits(b)
    api.lib.mm_b200_free_batch(b)
    one = api.opt_with(0)
    reads1, reads2 = _read_fq(r1), _read_fq(r2)
    assert len(got) == 2 * len(reads1)
    n_hits = 0
    for k in range(0, len(reads1), every):
        (n1, s1, _), (n2, s2, _) = reads1[k], reads2[k]
        want1, rep1 = api.map_frag(n1, [s1], one)
        want2, rep2 = api.map_frag(n2, [L.revcomp(s2) if flip2 else s2], one, len(s2) if flip2 else None)
        assert got[2 * k] == (want1[0], rep1), f"pair {k} mate 1"
        assert got[2 * k + 1] == (want2[0], rep2), f"pair {k} mate 2"
        n_hits += len(want1[0]) + len(want2[0])
    assert all(h[-1] == 0 for hits, _ in got for h in hits), "a hit has proper_frag set"
    return got, n_hits, list(pc)


@pytest.fixture(scope="module")
def synth(tmp_path_factory):
    if not (os.path.exists(SYN) and os.path.exists(NEW)):
        pytest.skip("needs build/mmsynth and build/minimap2-b200")
    d = tmp_path_factory.mktemp("nopair")
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "3000000", "3", "42"])
    subprocess.check_call([SYN, "sr", str(d / "ref.fa"), str(d / "r1.fq"), str(d / "r2.fq"), "4000", "46", "0.05"])
    _write_rc(d / "r2.fq", d / "r2rc.fq")
    return d


def test_api_sr_device_path(synth):
    api = Api(synth / "ref.fa", b"sr")
    try:
        got, n_hits, _ = _check_independent(api, synth / "r1.fq", synth / "r2.fq", True, every=4)
        assert n_hits > 1500
        # mm_b200_map_batches: several mini-batches, two in flight, each staged while the one before is mapped
        opt = api.opt_with(MM_F_INDEPEND_SEG)
        arr = (C.c_char_p * 2)(str(synth / "r1.fq").encode(), str(synth / "r2.fq").encode())
        reader = api.lib.mm_b200_open_reads(2, arr)
        bs = []
        while True:
            b = api.lib.mm_b200_read_batch(reader, C.byref(opt), 150_000)
            if not b:
                break
            bs.append(b)
        api.lib.mm_b200_close_reads(reader)
        assert len(bs) >= 6
        assert api.lib.mm_b200_map_batches(api.mi, C.byref(opt), 8, (C.c_void_p * len(bs))(*bs), len(bs), 0) == 0
        assert [x for b in bs for x in api.batch_hits(b)] == got
        for b in bs:
            api.lib.mm_b200_free_batch(b)
        # the joint mapping of the same pairs does pair them: the flag is what changed
        opt = api.opt_with(0)
        b = api.read_batch([synth / "r1.fq", synth / "r2.fq"], opt)
        assert api.lib.mm_b200_map_batch(api.mi, C.byref(opt), 8, b, 0) == 0
        joint = api.batch_hits(b)
        api.lib.mm_b200_free_batch(b)
        assert sum(h[-1] for hits, _ in joint for h in hits) > 1000
    finally:
        api.close()


def test_api_sr_paths_fixture(data):  # noqa: F811
    """re-chaining, warp hit trees, the heap replay and z-drop cuts under the flag: every pair is checked against the batch
    single-end path on r1 and revcomp(r2) (the same single-segment mapping as mm_map_frag, which checks every 8th pair)"""
    _write_rc(data / "r2.fq", data / "r2rc_np.fq")
    api = Api(data / "ref.fa", b"sr")
    try:
        L_ = api.lib
        got, n_hits, paths = _check_independent(api, data / "r1.fq", data / "r2.fq", True, every=8)
        assert n_hits > 1000
        one = api.opt_with(0)
        for fn, j in ((data / "r1.fq", 0), (data / "r2rc_np.fq", 1)):
            b = api.read_batch([fn], one)
            assert L_.mm_b200_map_batch(api.mi, C.byref(one), 8, b, 0) == 0
            want = api.batch_hits(b)
            L_.mm_b200_free_batch(b)
            reads = _read_fq(fn)
            for k, (w_hits, w_rep) in enumerate(want):
                if j == 1:  # back to the orientation of the read as it was read
                    ql = len(reads[k][1])
                    w_hits = [h[:3] + (ql - h[4], ql - h[3], 1 - h[5]) + h[6:] for h in w_hits]
                assert got[2 * k + j] == (w_hits, w_rep), f"pair {k} mate {j + 1}"
        # the batch under the flag: [0] rechained, [1] + [2] heap replays, [3] warp_tree, [4] zdrop_rounds, [5] zdrop_cuts.  Equal
        # positions in the seed merge come mostly from overlapping mates of one fragment, so the heap replay is rare here
        assert paths[0] > 100 and paths[3] > 100, paths
        assert paths[1] + paths[2] >= 1, paths
        assert paths[5] > 10 and paths[4] >= 1, paths
    finally:
        api.close()


def test_api_long_read_host_path(tmp_path):
    """-x map-ont --frag=yes on two files: the host stages (stage_hits / stage_finish); pe_ori = 0 flips nothing"""
    if not os.path.exists(SYN):
        pytest.skip("needs build/mmsynth")
    d = tmp_path
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "3000000", "3", "42"])
    subprocess.check_call([SYN, "long", str(d / "ref.fa"), str(d / "long.fq"), "120", "47", "4000"])
    reads = _read_fq(d / "long.fq")
    with open(d / "l1.fq", "wb") as f1, open(d / "l2.fq", "wb") as f2:
        for k in range(0, len(reads) - 1, 2):
            f1.write(_fastq(b"lp%d/1" % k, reads[k][1], reads[k][2]))
            f2.write(_fastq(b"lp%d/2" % k, reads[k + 1][1], reads[k + 1][2]))
    api = Api(d / "ref.fa", b"map-ont")
    try:
        api.opt.flag |= MM_F_FRAG_MODE
        assert api.opt.pe_ori == 0
        _, n_hits, _ = _check_independent(api, d / "l1.fq", d / "l2.fq", False)
        assert n_hits > 50
    finally:
        api.close()


def test_mm_map_frag_ignores_flag(synth):
    """the reference's mm_map_frag maps the segments it is given jointly whatever MM_F_INDEPEND_SEG says"""
    api = Api(synth / "ref.fa", b"sr")
    try:
        joint, indep = api.opt_with(0), api.opt_with(MM_F_INDEPEND_SEG)
        r1, r2 = _read_fq(synth / "r1.fq"), _read_fq(synth / "r2.fq")
        n_proper = 0
        for k in range(0, len(r1), 20):
            segs = [r1[k][1], L.revcomp(r2[k][1])]
            a = api.map_frag(r1[k][0], segs, joint)
            b = api.map_frag(r1[k][0], segs, indep)
            assert a == b, f"pair {k}"
            n_proper += sum(h[-1] for hits in a[0] for h in hits)
        assert n_proper > 50
    finally:
        api.close()


# ---------------------------------------------------------------------------------------------------- CLI

def _run(args, cwd):
    p = subprocess.run([NEW] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    return [l for l in p.stdout.decode().split("\n") if l and not l.startswith("@")]


def _by_read(lines):
    """records grouped by read, in order (each read's records are consecutive)"""
    out = []
    for l in lines:
        n = l.split("\t", 1)[0]
        if out and out[-1][0] == n:
            out[-1][1].append(l)
        else:
            out.append((n, [l]))
    return out


_PAIR_BITS = 0x1 | 0x2 | 0x8 | 0x20 | 0x40 | 0x80


def _toggle_sa(v):
    """SA:Z: value with every strand toggled"""
    out = []
    for e in v.split(";"):
        if e:
            x = e.split(",")
            x[2] = "+-"[x[2] == "+"]
            e = ",".join(x)
        out.append(e)
    return ";".join(out)


def _sam_norm(line, mate2):
    """a SAM record without its pairing fields; a mate-2 record of the paired run is brought to the single-end run on revcomp(r2)"""
    f = line.split("\t")
    name = f[0][:-2] if f[0][-2:] in ("/1", "/2") else f[0]
    flag = int(f[1]) & ~_PAIR_BITS
    if flag & 0x4:
        f[2], f[3] = "*", "0"  # an unmapped read is placed at its mate's primary in a pair
    if mate2:
        if not flag & 0x4:
            flag ^= 0x10
            for i in range(11, len(f)):
                if f[i].startswith("SA:Z:"):
                    f[i] = "SA:Z:" + _toggle_sa(f[i][5:])
        elif f[9] != "*":
            f[9] = L.revcomp(f[9].encode()).decode()
            f[10] = f[10][::-1]
    return "\t".join([name, str(flag)] + f[2:6] + f[9:])


def _paf_norm(line, l_seq=None):
    """a PAF record of the single-end run on revcomp(r2) in the read's own orientation (l_seq given), or as it is"""
    f = line.split("\t")
    if l_seq is not None:
        qs, qe = int(f[2]), int(f[3])
        f[2], f[3], f[4] = str(l_seq - qe), str(l_seq - qs), "+-"[f[4] == "+"]
    return "\t".join(f)


@pytest.mark.parametrize("extra", [[], ["--secondary=yes"], ["--cs", "--MD"], ["--paf"]], ids=lambda a: " ".join(a) or "sam")
def test_cli_equals_single_end(synth, extra):
    paf = extra == ["--paf"]
    x = ["-cx" if paf else "-ax", "sr"] + ([] if paf else extra) + ["-t", "8", "ref.fa"]
    got = _run(x[:2] + ["--no-pairing"] + x[2:] + ["r1.fq", "r2.fq"], synth)
    one1, one2 = _by_read(_run(x + ["r1.fq"], synth)), _by_read(_run(x + ["r2rc.fq"], synth))
    if paf:  # reads without a hit print nothing: pair the records by name
        d1, d2 = dict(one1), dict(one2)
        want = []
        for (n1, _, _), (n2, s2, _) in zip(_read_fq(synth / "r1.fq"), _read_fq(synth / "r2.fq")):
            want += d1.get(n1.decode(), []) + [_paf_norm(l, len(s2)) for l in d2.get(n2.decode(), [])]
        assert len(want) > 6000 and got == want
    else:
        assert len(one1) == len(one2) and len(one1) > 3000
        by = _by_read(got)  # paired QNAMEs are trimmed: a pair's records share one name
        assert len(by) == len(one1)
        for k, ((_, recs), (_, a), (_, b)) in enumerate(zip(by, one1, one2)):
            m1 = [_sam_norm(l, False) for l in recs if int(l.split("\t")[1]) & 0x40]
            m2 = [_sam_norm(l, True) for l in recs if int(l.split("\t")[1]) & 0x80]
            assert m1 == [_sam_norm(l, False) for l in a], f"pair {k} mate 1"
            assert m2 == [_sam_norm(l, False) for l in b], f"pair {k} mate 2"
            assert not any(int(l.split("\t")[1]) & 0x2 for l in recs)
    key = " ".join(["--no-pairing"] + x + ["r1.fq", "r2.fq"])
    if L.have_ref_bin():
        p = subprocess.run([L.REF_BIN_B] + x[:2] + ["--no-pairing"] + x[2:] + ["r1.fq", "r2.fq"], cwd=synth, stdout=subprocess.PIPE)
        assert p.returncode == 0
        want = [l for l in p.stdout.decode().split("\n") if l and not l.startswith("@")]
        assert len(want) == len(got)
        for i, (a, b) in enumerate(zip(want, got)):
            assert a == b, f"line {i}:\nref: {a[:300]}\nnew: {b[:300]}"
        return
    blob = "\n".join(got).encode()
    digest = {"bytes": len(blob), "sha256": hashlib.sha256(blob).hexdigest()}
    assert CLI_DIGESTS.get(key) == digest, f"{key!r}: {digest}"


def test_cli_two_gpus_same_bytes(synth):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    args = ["-ax", "sr", "--no-pairing", "-t", "8", "-K", "200k", "ref.fa", "r1.fq", "r2.fq"]
    assert _run(["--gpus", "2"] + args, synth) == _run(["--gpus", "1"] + args, synth)
