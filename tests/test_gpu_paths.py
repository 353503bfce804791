"""The kernels and code paths that only run for particular data must (a) actually run in the test suite and (b) give the
reference's bytes there.  The fixture is built for that: a 3 000-copy repeat family (minimizers between the two occurrence
cut-offs -> re-chain pass with thousands of chains per fragment), overlapping mates (equal positions meet in the seed merge),
reads with a block of mismatches (z-drop cuts), reads whose head is unrelated sequence (extension windows wider than the DP
band), and kilobase reads with an internal duplication mapped with the short-read preset (more merge lists than the rank
replay packs).  After each run the CLI's path counters / per-kernel launch counts (MM2_B200_PROFILE=1) are checked next to
the byte-for-byte comparison with oracle/_ref/minimap2_B, or with the output's digest recorded in tests/golden/digests.json where
the reference fork is not built."""
import os
import re
import subprocess
import numpy as np
import pytest
import _libs as L

pytestmark = pytest.mark.gpu
NEW = os.path.join(L.ROOT, "build", "minimap2-b200")


def _fastq(name, seq):
    return b"@" + name + b"\n" + seq + b"\n+\n" + b"I" * len(seq) + b"\n"


@pytest.fixture(scope="module")
def data(tmp_path_factory):
    if not os.path.exists(NEW):
        pytest.skip("needs build/minimap2-b200")
    d = tmp_path_factory.mktemp("paths")
    rng = np.random.default_rng(2024)
    ctg = [bytearray(L.rand_seq(rng, 2_000_000)) for _ in range(3)]
    elem = L.rand_seq(rng, 350)
    copies = []
    for i in range(3000):  # the high-copy family: every copy with its own 0-3 % divergence
        c, o = int(rng.integers(0, 3)), int(rng.integers(2000, 1_997_000))
        e = np.frombuffer(elem, dtype=np.uint8).copy()
        mut = rng.random(350) < rng.random() * 0.03
        e[mut] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, int(mut.sum()))]
        ctg[c][o:o + 350] = e.tobytes()
        copies.append((c, o))
    ctg = [bytes(c) for c in ctg]
    with open(d / "ref.fa", "wb") as f:
        for i, c in enumerate(ctg):
            f.write(b">chr%d\n" % (i + 1))
            f.write(b"\n".join(c[j:j + 80] for j in range(0, len(c), 80)) + b"\n")
    tr = bytes.maketrans(b"ACGT", b"CATG")
    r1, r2 = [], []

    def pair(name, frag, kind):
        if rng.random() < 0.5:
            frag = L.revcomp(frag)
        m1, m2 = bytearray(L.mutate(rng, frag[:150], 0.01, 0.0015, 0.0005)), bytearray(L.mutate(rng, L.revcomp(frag)[:150], 0.01, 0.0015, 0.0005))
        if kind == "zdrop" and len(m1) > 140:
            lo, ln = int(rng.integers(40, 70)), int(rng.integers(14, 45))
            m1[lo:lo + ln] = bytes(m1[lo:lo + ln]).translate(tr)
        if kind == "head" and len(m2) > 140:
            m2[:95] = L.rand_seq(rng, 95)
        r1.append(_fastq(name + b"/1", bytes(m1)))
        r2.append(_fastq(name + b"/2", bytes(m2)))

    for i in range(1200):  # fragments over a copy of the family
        c, o = copies[int(rng.integers(0, len(copies)))]
        st = o - int(rng.integers(20, 120))
        pair(b"rep%d" % i, ctg[c][st:st + int(rng.integers(300, 520))], "rep")
    for i in range(2500):  # unique sequence, short inserts: overlapping mates
        c = int(rng.integers(0, 3)); ins = int(np.clip(rng.normal(300, 70), 160, 600)); o = int(rng.integers(0, 2_000_000 - ins))
        pair(b"uni%d" % i, ctg[c][o:o + ins], ["uni", "uni", "uni", "zdrop", "head"][i % 5])
    open(d / "r1.fq", "wb").write(b"".join(r1))
    open(d / "r2.fq", "wb").write(b"".join(r2))
    with open(d / "kb.fq", "wb") as f:  # kilobase reads with an internal duplication, for the short-read preset single-end
        for i in range(24):
            c = int(rng.integers(0, 3)); o = int(rng.integers(0, 1_990_000))
            s = ctg[c][o:o + 2600]
            s = s[:1800] + s[600:1400] + s[1800:]
            f.write(_fastq(b"kb%d" % i, L.mutate(rng, s, 0.005, 0.001, 0.001)))
    with open(d / "long.fq", "wb") as f:
        for i in range(60):
            c = int(rng.integers(0, 3)); ln = int(rng.integers(1500, 9000)); o = int(rng.integers(0, 2_000_000 - ln))
            s = ctg[c][o:o + ln]
            f.write(_fastq(b"long%d" % i, L.mutate(rng, s if i % 2 else L.revcomp(s), 0.03, 0.03, 0.03)))
    return d


def _run(binary, args, cwd, profile=False):
    env = dict(os.environ, MM2_B200_PROFILE="1") if profile else None
    p = subprocess.run([binary] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    return [l for l in p.stdout.decode().split("\n") if not l.startswith("@PG")], p.stderr.decode()


def _stats(err):
    kern = {m.group(1): int(m.group(2)) for m in re.finditer(r"\[M::b200\] kernel (\S+)\s+(\d+) launches", err)}
    m = re.search(r"\[M::b200\] paths: (.*)", err)
    paths = {k: int(v) for k, v in re.findall(r"(\w+) (\d+)", m.group(1))} if m else {}
    return kern, paths


def _same_as_reference(args, got, cwd):
    if not L.have_ref_bin():
        L.check_digest("paths " + " ".join(args), got)
        return
    want, _ = _run(L.REF_BIN_B, args, cwd)
    assert len(want) == len(got)
    for i, (a, b) in enumerate(zip(want, got)):
        assert a == b, f"line {i}:\nref: {a[:300]}\nnew: {b[:300]}"
    L.record_reference_digest("paths " + " ".join(args), want)


def test_repeat_family_pairs(data):
    args = ["-ax", "sr", "-t", "8", "ref.fa", "r1.fq", "r2.fq"]
    got, err = _run(NEW, args, data, profile=True)
    _same_as_reference(args, got, data)
    kern, paths = _stats(err)
    assert paths.get("rechained", 0) > 100, paths            # the max_occ pass (map.c:353-375) and its CTA-per-fragment chain tail
    assert kern.get("k_chain_tail_block", 0) >= 1, kern
    assert paths.get("warp_tree", 0) > 100, paths             # hit trees of fragments with more than 32 chains
    assert paths.get("heap_rank_replay", 0) > 100, paths      # equal positions in the seed merge
    assert paths.get("zdrop_cuts", 0) > 10 and paths.get("zdrop_rounds", 0) >= 1, paths
    assert kern.get("k_ksw_tpj", 0) >= 1 and kern.get("k_ksw_dpx", 0) >= 1, kern   # both DP forms


def test_kilobase_reads_short_read_preset(data):
    args = ["-ax", "sr", "-t", "4", "ref.fa", "kb.fq"]
    got, err = _run(NEW, args, data, profile=True)
    _same_as_reference(args, got, data)
    kern, paths = _stats(err)
    assert paths.get("heap_literal_replay", 0) + paths.get("heap_rank_replay", 0) >= 1, paths


def test_long_reads_wavefront_dp(data):
    args = ["-ax", "map-ont", "-t", "8", "ref.fa", "long.fq"]
    got, err = _run(NEW, args, data, profile=True)
    _same_as_reference(args, got, data)
    kern, _ = _stats(err)
    assert kern.get("k_ksw_wave", 0) >= 1, kern
